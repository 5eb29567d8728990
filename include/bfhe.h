/*
 * bfhe.h -- C ABI of the B200-native gate-bootstrapping engine.
 *
 * This is the drop-in boundary beneath the reference's circuit evaluator.  Each entry point
 * names the lbcrypto::BinFHEContext call (and the call site in /root/reference) it replaces.
 * Plain pointers and sizes only; no C++ or torch types.  All functions return 0 on success and
 * a negative code on error (text from bfhe_last_error()); nothing throws across this boundary.
 *
 * Ciphertexts: an LWE ciphertext mod q is ct_words = n+1 uint32 words (a_0..a_{n-1}, b) stored in a
 * row of ct_stride words (ct_words rounded up to a multiple of 4).  A "slab" is a device array of
 * such rows; gates name their operands by row index, exactly like the reference's registers
 * (R<k> in the .out format, src/circuit.cpp:144-294).
 *
 * There is NO CPU fallback: every Eval* entry point runs hand-written sm_100a kernels and fails
 * with BFHE_ERR_CUDA when no device is available.
 */
#ifndef BFHE_H
#define BFHE_H
#include <stddef.h>
#include <stdint.h>
#ifdef __cplusplus
extern "C" {
#endif

/* enum values follow OpenFHE 1.0.x binfhe-constants.h (lbcrypto::BINFHE_PARAMSET / BINFHE_METHOD / BINGATE);
 * the reference only ever passes TOY / STD128_OPT and AP / GINX (src/circuit.cpp:69-86, src/utils.cpp:165-190) */
enum { BFHE_TOY = 0, BFHE_STD128_OPT = 5 };
enum { BFHE_AP = 0, BFHE_GINX = 1 };
enum { BFHE_OR = 0, BFHE_AND = 1, BFHE_NOR = 2, BFHE_NAND = 3, BFHE_XOR_FAST = 4, BFHE_XNOR_FAST = 5,
       BFHE_XOR = 6, BFHE_XNOR = 7, /* composite OR(AND(a,!b),AND(!a,b)) as src/gate.cpp:198-202 */
       BFHE_BOOTSTRAP = 8 /* BinFHEContext::Bootstrap: in1 ignored */ };
#define BFHE_NEG0 0x100u /* operand 0 passes through EvalNOT first (fused, no bootstrap) */
#define BFHE_NEG1 0x200u

enum { BFHE_OK = 0, BFHE_ERR_ARG = -1, BFHE_ERR_STATE = -2, BFHE_ERR_CUDA = -3, BFHE_ERR_FORMAT = -4,
       BFHE_ERR_ALIAS = -5 /* EvalBinGate(ct, ct): OpenFHE throws, src/gate.cpp:134 catches */,
       BFHE_ERR_NCCL = -6, BFHE_ERR_IO = -7 };

typedef struct {
  uint32_t paramset, method;
  uint32_t n, N, q;
  uint64_t Q, qKS;
  uint32_t baseKS, dKS, baseG, dG, baseR, dR;
  uint32_t ct_words, ct_stride;
} bfhe_params;

/* one gate of a wavefront: replaces one Gate::Evaluate task (src/gate.cpp:49, src/circuit.cpp:698-710) */
typedef struct {
  uint32_t op; /* BFHE_<gate> | BFHE_NEG0 | BFHE_NEG1 */
  uint32_t in0, in1, out; /* slab rows */
} bfhe_gate;

typedef struct bfhe_ctx bfhe_ctx;

/* ---- context: BinFHEContext::GenerateBinFHEContext(set, method)  (src/circuit.cpp:88) ---- */
bfhe_ctx *bfhe_create(int paramset, int method, int device /* CUDA ordinal, -1 = host-only (keygen/encrypt/decrypt) */);
void bfhe_destroy(bfhe_ctx *);
int bfhe_get_params(const bfhe_ctx *, bfhe_params *out);
const char *bfhe_last_error(void);
/* launch stream for every subsequent kernel: a cudaStream_t (e.g. torch's current stream; NULL = the legacy default
 * stream), or use_own != 0 to go back to the context's private non-blocking stream (the initial state) */
int bfhe_set_stream(bfhe_ctx *, void *cuda_stream, int use_own);
int bfhe_sync(bfhe_ctx *);

/* ---- keys: KeyGen() / BTKeyGen(sk)  (src/circuit.cpp:90-91) ----
 * Randomness contract (keygen, btkeygen, encrypt, circuit_set_input): every secret, mask and noise term is drawn from a ChaCha20
 * stream.  seed == 0 keys the stream with 256 bits of OS entropy (getrandom): the secure default, equivalent to OpenFHE's self-seeding
 * PRNG that the reference relies on.  seed != 0 derives the stream from the 64-bit seed alone: reproducible keys / ciphertexts for
 * tests, oracle parity and benchmarks, and therefore NOT confidential.  For sharded (multi-rank) evaluation generate the keys on one
 * rank with seed 0 and distribute the blob (bfhe_export_keys -> broadcast -> bfhe_import_keys); do not share a constant seed. */
int bfhe_keygen(bfhe_ctx *, uint64_t seed);   /* LWE secret key (host) */
int bfhe_btkeygen(bfhe_ctx *, uint64_t seed); /* bootstrapping + key-switching keys (host), uploaded if a device is attached */
/* flat key blob ("same serialized keys" contract, SURVEY 5 checkpoint/resume): layout documented in DESIGN.md:
 *   header{magic "BFHEKEY1", version, params, has_sk, ksk_elem_bytes, Q, qKS, bk_words, ksk_elems}
 *   sk[n] int32 | BK coefficient form uint32 | KSK [N][baseKS][dKS][n+1] uint16 (qKS<=2^16) or uint32 */
size_t bfhe_keyblob_size(const bfhe_ctx *);
int bfhe_export_keys(const bfhe_ctx *, void *buf, size_t cap, int include_sk);
/* either blob, BFHEKEY1 or BFHEKEY2 (below); the parameters must match this context, else BFHE_ERR_FORMAT */
int bfhe_import_keys(bfhe_ctx *, const void *buf, size_t len);
int bfhe_save_keys(const bfhe_ctx *, const char *path, int include_sk);
int bfhe_load_keys(bfhe_ctx *, const char *path);

/* ---- compact evaluation keys: the public masks come from a seed ----
 * Most of a key blob is uniform masks that carry no secret: n of the n+1 words of every KSK row, and column 0 of every RGSW row of the
 * BK.  bfhe_btkeygen_compact generates the same kinds of keys as bfhe_btkeygen, with the same noise, and leaves the context in the same
 * state, but every mask is the expansion of a 256-bit public MASK SEED that the context keeps.  Its blob, BFHEKEY2, then carries only the
 * seed and the bodies: at STD128_OPT about 33.4 MB instead of 329.5 MB (GINX) and 1.02 GB instead of 2.30 GB (AP).
 *   mask seed: seed == 0 -> 256 bits of OS entropy, drawn independently of the secret stream; seed != 0 -> 256 bits of a dedicated stream
 *              of the secret SeedKey (reproducible for tests, and ChaCha20 output reveals nothing about its key).
 *   expansion: mask row r is the ChaCha20 keystream (RFC 8439 block function, 64-bit block counter from 0 in words 12-13, 64-bit nonce
 *              in words 14-15) with key = mask seed (eight little-endian words) and nonce = r.  Coefficient t of the row is the
 *              little-endian 128-bit integer of keystream words 4t .. 4t+3, reduced mod the row's modulus m (qKS for the KSK, Q for the
 *              BK): statistical distance from uniform below m / 2^128 per coefficient, no rejection, so one ChaCha block gives four
 *              coefficients and any of them can be computed alone.
 *   rows:      KSK row (i, j, k) (i < N, digit value j < baseKS, digit k < dKS) is r = (i * baseKS + j) * dKS + k; BK mask polynomial p is
 *              r = 2^40 + p, where p counts the column-0 polynomials in BFHEKEY1 order (RGSW t, row l: p = t * 2dG + l).
 *   bodies:    KSK b = <a,s> + e + z_i * j * baseKS^k mod qKS, as bfhe_btkeygen.  BK row l of an RGSW of m (m = 1 or 0 for GINX,
 *              +-X^mm for AP): odd rows b = a*z + e + m*g^(l/2), as bfhe_btkeygen; even rows, whose message bfhe_btkeygen adds to the
 *              mask, b = a*z + e - m*g^(l/2)*z, so the public mask never carries the message.  The phase b - a*z is unchanged, and the
 *              kernels see an ordinary RGSW key.
 * SECURITY: the mask seed is public.  It is drawn fresh by every call, so two key sets never share one; never reuse a mask seed for
 * another key set (two key sets with one seed and different secrets would share their masks).
 * Layout of BFHEKEY2: the BFHEKEY1 header with magic "BFHEKEY2", version 1 (the same fields and values) | mask seed, 32 bytes |
 *   sk[n] int32 (zero without the secret key) | BK bodies: the column-1 polynomials in BFHEKEY1 order, coefficient form, uint32 |
 *   KSK bodies [N][baseKS][dKS], uint16 when qKS <= 2^16 else uint32; each section padded to 8 bytes, as in BFHEKEY1.
 * Import checks every body word against its modulus (BFHE_ERR_FORMAT naming the section and index, before any device work, leaving the
 * previous keys in place).  A device context uploads the bodies and generates the masks on the GPU; it keeps the bodies, not the full
 * keys, on the host, and bfhe_export_keys / bfhe_export_openfhe_json expand them on the host when called.  A host-only context expands
 * them on import. */
int bfhe_btkeygen_compact(bfhe_ctx *, uint64_t seed);
size_t bfhe_keyblob_compact_size(const bfhe_ctx *);
/* BFHE_ERR_STATE when the keys have no mask seed (bfhe_btkeygen, a BFHEKEY1 import, an OpenFHE JSON import) */
int bfhe_export_keys_compact(const bfhe_ctx *, void *buf, size_t cap, int include_sk);

/* ---- compact fresh ciphertexts: a client's inputs as a public mask seed and one body word per bit ----
 * n of the n+1 words of a fresh encryption are its uniform mask, which carries no secret.  bfhe_encrypt_compact draws every mask from a
 * public seed, so the blob, BFHECTS1, holds that seed and one body per bit: an AES-128 block (256 bits) is 576 bytes instead of 516 KB of
 * full rows at STD128_OPT.  Only fresh encryptions can be compact; bootstrapped ciphertexts and the evaluator's outputs stay full rows.
 *   mask seed: 256 bits, fresh on every call.  seed == 0 -> OS entropy, independent of the secret stream; seed != 0 -> a dedicated stream
 *              of the secret SeedKey (reproducible and not confidential, as for every nonzero seed; a different stream from the mask
 *              seed of bfhe_btkeygen_compact).
 *   expansion: row g (g = 0 .. count-1) has mask row r = g under this seed, by the rule of the compact keys above: ChaCha20 keyed with the
 *              seed, nonce r, coefficient t = keystream words 4t .. 4t+3 as a little-endian 128-bit integer mod q.  q is a power of two,
 *              so the reduction is exact and uniform.
 *   body:      b_g = <a_g, s> + e_g + (bits[g] % 4) * q/4 mod q, the message convention of bfhe_encrypt; e_g is the Gaussian noise of
 *              bfhe_encrypt drawn from stream 2^48 + g of the secret SeedKey (a range no other call uses).
 * Layout of BFHECTS1, little-endian: 64-byte header {magic "BFHECTS1", u32 version = 1, u32 paramset, u32 n, u32 q, u64 count, the 32-byte
 *   mask seed} | count uint16 bodies, zero-padded to 8 bytes.  Size 64 + pad8(2 * count).
 * Every reader checks on the host, before any device work, and answers BFHE_ERR_FORMAT naming what failed: magic and version; paramset,
 *   n and q equal to the context's; the exact length; every body below q (naming the first bad index); zero padding bytes.
 * SECURITY: the mask seed is public and the noise comes only from the secret stream.  Never reuse a mask seed for a second batch under
 * the same key: identical masks expose the differences of the messages.  bfhe_encrypt_compact draws a new one on every call. */
size_t bfhe_ct_compact_size(const bfhe_ctx *, size_t count);
/* on the host, with the secret key (BFHE_ERR_STATE without it); works on host-only contexts.  blob holds bfhe_ct_compact_size bytes. */
int bfhe_encrypt_compact(const bfhe_ctx *, const uint8_t *bits, size_t count, uint64_t seed, void *blob, size_t cap);
/* the blob's count full rows of ct_stride words (padding words zero) into cts (cap_rows rows).  on_device == 0: host memory, works on any
 * context, with or without keys.  on_device != 0: memory of the context's device, 16-byte aligned (else BFHE_ERR_ARG), written by one
 * expansion launch on the launch stream; returns after the rows are written.  A host-only context gives BFHE_ERR_CUDA. */
int bfhe_expand_cts(bfhe_ctx *, const void *blob, size_t len, uint32_t *cts, size_t cap_rows, int on_device);

/* ---- OpenFHE 1.0.x object exchange (SURVEY 8 row f-3; the reference's crypto is find_package(OpenFHE), CMakeLists.txt:8, "Tested with
 * OpenFHE v.1.0.1", Release_Notes.md:4) ----
 * cereal JSON archives as OpenFHE's own Serial::SerializeToFile(path, obj, SerType::JSON) writes them (the reference itself never
 * serialises): the LWE secret key (LWEPrivateKey), the refresh key (cc.GetRefreshKey(), RingGSWACCKey), the switching key
 * (cc.GetSwitchKey(), LWESwitchingKey) and single LWE ciphertexts.  Refresh-key polynomials are taken in EVALUATION format (OpenFHE's
 * order: Cooley-Tukey bit-reversed, smallest primitive 2N-th root) or COEFFICIENT format, per polynomial as its "f" member says.
 * Importing both the refresh and the switching key leaves the context exactly as after bfhe_btkeygen.  A file whose ring modulus is
 * not this context's Q is refused with BFHE_ERR_FORMAT (DESIGN.md section 3).  The layout is restated from the 1.0.x sources from
 * memory -- OpenFHE is not available in this build environment -- so parity against a real OpenFHE file is UNPINNED until a
 * maintainer runs tools/openfhe_export_keys.cpp (INTEGRATION.md "Closing the parity gap").  cereal's portable-binary form is
 * positional and cannot be checked offline; it is deliberately not offered. */
enum { BFHE_OFHE_SECRET_KEY = 0, BFHE_OFHE_REFRESH_KEY = 1, BFHE_OFHE_SWITCH_KEY = 2 };
int bfhe_import_openfhe_json(bfhe_ctx *, int what, const char *path);
int bfhe_export_openfhe_json(const bfhe_ctx *, int what, const char *path);
int bfhe_import_openfhe_ct_json(const bfhe_ctx *, const char *path, uint32_t *ct_row /* ct_stride words */);
int bfhe_export_openfhe_ct_json(const bfhe_ctx *, const uint32_t *ct_row, const char *path);

/* ---- host-side LWE: Encrypt(sk, bit, FRESH) / Decrypt(sk, ct, &res)  (src/circuit.cpp:506,800; src/gate.cpp:72..) ---- */
int bfhe_encrypt(const bfhe_ctx *, const uint8_t *bits, size_t count, uint64_t seed, uint32_t *ct_host /* count*ct_stride */);
int bfhe_decrypt(const bfhe_ctx *, const uint32_t *ct_host, size_t count, uint8_t *out /* floor(4r/q) in 0..3 */);

/* ---- device slabs (wire storage; replaces Wire::ct shared_ptrs, src/wire.h:46-73) ---- */
int bfhe_slab_alloc(bfhe_ctx *, size_t rows, uint32_t **dev_ptr);
int bfhe_slab_free(bfhe_ctx *, uint32_t *dev_ptr);
int bfhe_slab_upload(bfhe_ctx *, uint32_t *dev_slab, size_t first_row, const uint32_t *host, size_t rows);
int bfhe_slab_download(bfhe_ctx *, const uint32_t *dev_slab, size_t first_row, uint32_t *host, size_t rows);

/* ---- the hot path ---- */
/* EvalNOT(ct) for a batch (src/gate.cpp:112) */
int bfhe_eval_not_batch(bfhe_ctx *, uint32_t *dev_slab, const uint32_t *in_rows, const uint32_t *out_rows, size_t count);
/* EvalBinGate(gate, ct1, ct2) for one wavefront of independent gates (src/gate.cpp:133,146,172,200-202).
 * gates is a HOST array; XOR/XNOR expand to the reference's 3-bootstrap composite.  Asynchronous on the stream. */
int bfhe_eval_bingate_batch(bfhe_ctx *, uint32_t *dev_slab, const bfhe_gate *gates, size_t count);
/* Bootstrap(ct) for a batch (what Encrypt's BOOTSTRAPPED default applies to every input, src/circuit.cpp:506) */
int bfhe_bootstrap_batch(bfhe_ctx *, uint32_t *dev_slab, const uint32_t *in_rows, const uint32_t *out_rows, size_t count);
/* end-to-end form with HOST buffers: H2D of the input slab rows, the wavefront, D2H of the produced rows.
 * in_host holds rows [0, in_rows) of the slab; gate.out rows are >= in_rows and < in_rows + out_rows.  The padding words of every
 * output row are zero.
 * Concurrent calls on one context may be combined into one wave: a call that finds no batch in flight launches at once with whatever
 * is queued; calls that arrive while a batch runs queue up and go together as the next batch.  Results are identical to separate calls
 * (a gate's words do not depend on the batch it ran in), and each call returns after its own rows are written.  Each call's arguments
 * (pointers, row ranges, op, the alias rule) are checked in its own thread before it joins, so a bad call fails alone; a CUDA failure
 * during a batch fails every call in it, each with the message in its own bfhe_last_error(). */
int bfhe_eval_bingate_host(bfhe_ctx *, const bfhe_gate *gates, size_t count, const uint32_t *in_host, size_t in_rows,
                           uint32_t *out_host, size_t out_rows);
/* EvalNOT(ct) on the host, for count rows of HOST memory: needs no device and works on host-only contexts.  The words of the device
 * EvalNOT: a_i -> (q - a_i) mod q, b -> (q/4 + q - b) mod q; padding words are written as zero.  Every input word a_0 .. a_{n-1}, b
 * must be below q, else BFHE_ERR_FORMAT naming the first bad row, and nothing is written.  ct_out may equal ct_in. */
int bfhe_eval_not_host(const bfhe_ctx *, const uint32_t *ct_in, size_t count, uint32_t *ct_out);

/* ---- measurement hooks ---- */
/* when enabled, every hot-path launch is bracketed by CUDA events on the launch stream */
int bfhe_profile_enable(bfhe_ctx *, int on);
/* kernel: 0 = blind rotation, 1 = key switch, 2 = EvalNOT; returns accumulated device ms and launch count, then resets */
int bfhe_profile_read(bfhe_ctx *, int kernel, double *ms, uint64_t *launches);
/* integer-pipe microbenchmark: measured 32-bit multiply-class instructions/s (IMAD, IMAD.HI, IMAD.WIDE) */
int bfhe_microbench_int(bfhe_ctx *, int which, double *ginstr_per_s);

/* ---- stage-level entry points (parity tests against the oracle; same kernels the hot path launches) ---- */
int bfhe_dbg_ntt_roundtrip(bfhe_ctx *, const uint32_t *poly_host, size_t npoly, uint32_t *fwd_inv_host, uint32_t *prod_host,
                           const uint32_t *poly2_host);
/* blind rotation only: acc in coefficient form (2N words per gate) */
int bfhe_dbg_blind_rotate(bfhe_ctx *, uint32_t *dev_slab, const bfhe_gate *gates, size_t count, uint32_t *acc_host);
/* test hook: force the blind-rotation form.  0 = cost model; 1, 2, 4 = that many gates per CTA (first-generation throughput
 * kernel); 8 = one gate per CTA, TMA-staged key (latency kernel); 32 = one gate on a 2-CTA thread-block cluster (STD128_OPT GINX);
 * 128 = one gate on a slot-sliced 4-CTA cluster (STD128_OPT, GINX and AP).  16 and 64 named round-1 forms that no longer exist. */
int bfhe_dbg_set_gates_per_cta(bfhe_ctx *, int gates_per_cta);
/* how many gates the 2-CTA / 4-CTA cluster forms keep co-resident on this device (cudaOccupancyMaxActiveClusters; differs between GPUs) */
int bfhe_dbg_cluster_limits(bfhe_ctx *, int *cl2_gates, int *cl4_gates);
/* imports a BFHEKEY2 blob as bfhe_import_keys does on a device context (same kernels and buffers) and writes the BFHEKEY1 blob the device
 * expansion produced: the BK staging buffer as downloaded, the device KSK restored to [N][baseKS][dKS][n+1] on the host.  full_blob holds
 * bfhe_keyblob_size bytes; the context keeps the imported keys. */
int bfhe_dbg_expand_keys(bfhe_ctx *, const void *compact_blob, size_t len, void *full_blob, size_t cap);
/* test hook for the combining of bfhe_eval_bingate_host: while hold != 0, calls queue and nothing launches, not even from an idle
 * context; hold = 0 launches everything queued as one batch (in one of the waiting callers' threads).  Returns the number of calls
 * that were queued when it was called (>= 0), so a test can wait until every caller has joined, or BFHE_ERR_ARG. */
int bfhe_dbg_hold_batches(bfhe_ctx *, int hold);

/* ---- circuit evaluator: mirrors class Circuit (src/circuit.h:56-72), level-synchronous ---- */
typedef struct bfhe_circuit bfhe_circuit;
bfhe_circuit *bfhe_circuit_create(bfhe_ctx *);
void bfhe_circuit_destroy(bfhe_circuit *);
int bfhe_circuit_read_file(bfhe_circuit *, const char *path);             /* Circuit::ReadFile (.out assembler format) */
int bfhe_circuit_read_bristol(bfhe_circuit *, const char *path, int new_format); /* analyze+assemble without the text round trip */
/* netlist from arrays / back to arrays / emitted as the reference's ".out" text.  kind[] uses GateEnum order
 * {INPUT, OUTPUT, NOT, AND, OR, XOR, DFF, LUT3, LUT4} (src/gate.h:51), then the native single-bootstrap gate types of EvalBinGate and
 * the composite XNOR: {NAND, NOR, XNOR, XOR_FAST, XNOR_FAST}.  INPUT: in0 = bus, in1 = bit, out = wire; OUTPUT: in0 = wire, out = bit;
 * DFF: in0 = D, out = Q (state 0 after Reset; Clock() may be called repeatedly, each call latches D -- the reason the reference's
 * method is called Clock(), README.md:55); LUT3 / LUT4 (stubs in the reference, src/gate.cpp:220-225): in0..in3 and a truth table whose
 * bit (in0 | in1 << 1 | in2 << 2 | in3 << 3) is the output, lowered at load to <= 5 / <= 13 two-input gates (_ex entry point).
 * ".out" grammar of the additions: "R3 = NAND(R1, R2)", "R5 = DFF(R4)", "R9 = LUT3(R1, R2, R3, 0xE8)", "R9 = LUT4(R1, R2, R3, R4, 0x6996)". */
int bfhe_circuit_load_netlist(bfhe_circuit *, const uint8_t *kind, const uint32_t *in0, const uint32_t *in1, const uint32_t *out,
                              size_t count, uint32_t n_wires, const uint32_t *in_bits, uint32_t n_in_buses, uint32_t out_bits);
int bfhe_circuit_load_netlist_ex(bfhe_circuit *, const uint8_t *kind, const uint32_t *in0, const uint32_t *in1, const uint32_t *in2,
                                 const uint32_t *in3, const uint32_t *table, const uint32_t *out, size_t count, uint32_t n_wires,
                                 const uint32_t *in_bits, uint32_t n_in_buses, uint32_t out_bits);
int bfhe_circuit_get_netlist(const bfhe_circuit *, uint8_t *kind, uint32_t *in0, uint32_t *in1, uint32_t *out, size_t cap,
                             uint32_t *count, uint32_t *n_wires);
int bfhe_circuit_write_out(const bfhe_circuit *, const char *path);
int bfhe_circuit_set_flags(bfhe_circuit *, int plaintext, int encrypted, int verify); /* setPlaintext/Encrypted/Verify */
int bfhe_circuit_info(const bfhe_circuit *, uint32_t *n_inputs, uint32_t *input_bits /*[8]*/, uint32_t *n_output_bits,
                      uint32_t *n_gates, uint32_t *n_bootstraps, uint32_t *n_levels, uint32_t *max_width);
/* multi-GPU: shard every level over world ranks; comm_id = 128-byte ncclUniqueId distributed by the caller.  From here on set_sharding,
 * set_wave_capacity, set_shard_threshold, set_flags, set_input and clock are COLLECTIVE: every rank makes the same calls in the same order
 * (they exchange launch costs and memory handles, and a rank's Clock stores into its peers' slabs) */
int bfhe_circuit_set_sharding(bfhe_circuit *, int rank, int world, const void *nccl_unique_id);
int bfhe_get_nccl_unique_id(void *out128);
/* how the ranks exchange a sharded level's output ciphertexts: 0 = single rank; 2 = the key-switch kernel stores every output into every
 * rank's slab itself (peer slabs mapped with CUDA IPC, stores over NVLink, one flag per rank and level -- chosen when every rank could
 * map every slab); 1 = one ncclAllGather per level (fallback, or BFHE_EXCHANGE=nccl in the environment).  Valid after the first
 * encrypted SetInput. */
int bfhe_circuit_exchange_mode(const bfhe_circuit *);
/* schedule: 0 = the reference's ASAP waves (src/circuit.cpp:593-677), one launch per level; n > 0 = ready gates packed into
 * waves of at most n bootstraps by longest remaining path; -1 (default) = one gate per SM and rank when a device is attached,
 * ASAP otherwise.  Ciphertexts do not depend on the schedule.  bfhe_circuit_info always reports the ASAP statistics. */
int bfhe_circuit_set_wave_capacity(bfhe_circuit *, int max_bootstraps_per_wave);
/* multi-GPU: levels with fewer than min_bootstraps bootstraps are computed redundantly by every rank and skip the exchange
 * (SURVEY 8(e)); 0 = shard every level; -1 (default) = per level by the measured cost model (device attached), else shard all */
int bfhe_circuit_set_shard_threshold(bfhe_circuit *, int min_bootstraps);
int bfhe_circuit_reset(bfhe_circuit *);                                     /* Circuit::Reset */
int bfhe_circuit_set_input(bfhe_circuit *, const uint8_t *bits, size_t nbits, uint64_t seed); /* Circuit::SetInput (all input buses concatenated) */
int bfhe_circuit_clock(bfhe_circuit *, uint8_t *out_bits, size_t cap, uint8_t *plain_out_bits); /* Circuit::Clock */
/* ---- evaluation with the evaluation keys only (a context that imported bfhe_export_keys(..., include_sk = 0)) ----
 * Circuit::SetInput on ciphertexts.  Needs evaluation keys only, never the secret key.  cts: nbits rows of ct_stride words, the input
 * buses concatenated in SetInput's bit order; on_device != 0: memory on the context's device, read in order on the launch stream
 * (bfhe_set_stream), else host memory.  Level 0 bootstraps them, exactly as it bootstraps SetInput's fresh encryptions.
 * Input contract: every word a_0 .. a_{n-1}, b is below q, else BFHE_ERR_FORMAT naming the first bad row, and the circuit is left
 * without input (Clock fails with BFHE_ERR_STATE until the next SetInput).  Padding words are ignored and stored as zero.
 * Modes: encrypted mode with plaintext and verify mode off, else BFHE_ERR_STATE (ciphertext inputs have no plaintext).  Argument and
 * state errors are reported before the device is touched.
 * Flip-flops power up from the trivial encryption of 0 (all-zero row), bootstrapped into the latch row: they decrypt exactly as after
 * SetInput(bits), whose power-up value is Encrypt(0), but the state rows' ciphertexts differ.
 * Sharded circuits (world > 1): collective; rank 0's rows are used and broadcast with rank 0's validation status, so every rank returns
 * the same code.  Other ranks may pass NULL.
 * After this call bfhe_circuit_clock (bits) decrypts as usual when the context holds the secret key, and fails with BFHE_ERR_STATE
 * before launching anything when it does not. */
int bfhe_circuit_set_input_ct(bfhe_circuit *, const uint32_t *cts, size_t nbits, int on_device);
/* bfhe_circuit_set_input_ct from a BFHECTS1 blob (bfhe_encrypt_compact): the masks are generated on the GPU straight into the circuit's
 * fresh input rows.  Modes, flip-flop power-up and the "without input on error" rule are those of bfhe_circuit_set_input_ct.  The blob's
 * checks give BFHE_ERR_FORMAT; count != the circuit's input bits gives BFHE_ERR_ARG.  Sharded circuits: collective; only rank 0's blob is
 * read (other ranks may pass NULL), and a blob rank 0 refuses still goes through the broadcast, so every rank returns the same code. */
int bfhe_circuit_set_input_compact(bfhe_circuit *, const void *blob, size_t len);
/* Circuit::Clock with the outputs left encrypted: out_bits rows of ct_stride words (padding words zero) into out_cts, host or device
 * memory (on_device as above).  An output that reads its wire through NOT comes out as EvalNOT of that row, so it decrypts to what
 * bfhe_circuit_clock returns.  Encrypted mode without verify mode; works after either SetInput form and needs no secret key.  Every rank
 * of a sharded circuit returns all outputs.  Returns after the rows are written. */
int bfhe_circuit_clock_ct(bfhe_circuit *, uint32_t *out_cts, size_t cap_rows, int on_device);
int bfhe_circuit_stats(const bfhe_circuit *, double *device_ms, double *host_ms, uint64_t *verify_mismatches);
/* the schedule in use: wave capacity (0 = ASAP), levels incl. the input-bootstrap level, levels that are sharded, and the four launch
 * costs (ms: 4-CTA cluster, 2-CTA cluster, one gate per SM, four gates per SM) the planner used -- measured by a start-up probe on the
 * first encrypted SetInput when the capacity is left to the cost model */
int bfhe_circuit_get_schedule(const bfhe_circuit *, uint32_t *wave_cap, uint32_t *n_levels, uint32_t *n_sharded, double *cost_ms4);
/* per-level plan, for tests of the sharding logic: gates of level L assigned to `rank` of `world`; *rows_per_rank == 0 with
 * world > 1 means the level is not sharded (every rank evaluates all of it, no exchange follows) */
int bfhe_circuit_level_plan(const bfhe_circuit *, uint32_t level, int rank, int world, bfhe_gate *out, size_t cap,
                            uint32_t *count, uint32_t *first_row, uint32_t *rows_per_rank);
/* plan internals for tests: total slab rows, first fresh-encryption row, level count incl. the input-bootstrap
 * level 0, slab row of every output bit (bit 31 set = read through NOT), and the EvalNOT pairs of one level */
int bfhe_circuit_plan_misc(const bfhe_circuit *, uint32_t *total_rows, uint32_t *fresh_base, uint32_t *n_levels_incl_input,
                           uint32_t *out_rows, uint32_t *not_count, uint32_t level, uint32_t *not_pairs);
int bfhe_circuit_use_graph(bfhe_circuit *, int on); /* one CUDA graph per circuit instead of per-level launches (default on) */
int bfhe_circuit_download_slab(bfhe_circuit *, uint32_t *host, size_t rows_cap); /* every wire ciphertext, for parity tests */
int bfhe_circuit_dump_gate_count(const bfhe_circuit *, uint32_t *in, uint32_t *out, uint32_t *and_, uint32_t *or_,
                                 uint32_t *xor_, uint32_t *not_);
int bfhe_circuit_dump_gate_count_ex(const bfhe_circuit *, uint32_t *counts8 /* DFF, LUT3, LUT4, NAND, NOR, XNOR, XOR_FAST, XNOR_FAST */);
/* Circuit::dumpNetList (what = 0: wire name -> names of the gates reading it, in the reference's map order) / Circuit::dumpGates
 * (what = 1: input gate names, then all gate names) as text (src/circuit.cpp:844-865); *needed = length without the final 0 */
int bfhe_circuit_dump_text(const bfhe_circuit *, int what, char *buf, size_t cap, size_t *needed);
/* clocked circuits, for tests of the plan: per flip-flop {row D is read from | bit 31 = through EvalNOT, state row (Q), latch row,
 * row of the fresh Encrypt(0) that the first clock after Reset bootstraps into the latch row} */
int bfhe_circuit_dff_plan(const bfhe_circuit *, uint32_t *n_dff, uint32_t *quads, size_t cap_dffs);

#ifdef __cplusplus
}
#endif
#endif
