--[[ ganrev.lua -- LuaJIT-FFI binding of libganrev_cuda.so (include/ganrev.h).

Drop-in arithmetic for aleju/gan-reverser's apply_r.lua: the models.lua G/R constructors and
apply_r.lua's search, cluster, fix and anomaly modes keep their names and call this module
instead of nn / cudnn / unsup / torch.dist.  No cutorch, no cudnn, no CPU fallback.

NOT EXECUTED IN THIS REPOSITORY'S CI: the build image has no lua/luajit/th.  Every call below
is mirrored one-to-one by gan-reverser_b200/_lib.py (ctypes), which is what the tests drive.

Usage (see INTEGRATION.md):
    local ganrev = require 'ganrev'
    local ctx = ganrev.new(OPT.gpu)                       -- replaces cutorch.setDevice(OPT.gpu + 1)
    MODEL_G = ganrev.wrap_G(ctx, tmp.G, {1, 32, 32}, 100)  -- flattens the trained nn.Sequential
    images  = MODEL_G:forward(noise)
]]
local ffi = require 'ffi'
require 'torch'

ffi.cdef[[
int usleep(unsigned int usec);
typedef struct ganrev_ctx ganrev_ctx;
int         ganrev_version(void);
int         ganrev_create(ganrev_ctx** out, int device);
void        ganrev_destroy(ganrev_ctx* ctx);
const char* ganrev_last_error(const ganrev_ctx* ctx);
int ganrev_comm_unique_id(ganrev_ctx* ctx, void* out, size_t cap, size_t* len);
int ganrev_comm_init(ganrev_ctx* ctx, int world, int rank, const void* uid, size_t len);
int ganrev_load_G(ganrev_ctx* ctx, int C, int H, int W, int noise_dim, const float* blob, size_t n_floats);
int ganrev_load_R(ganrev_ctx* ctx, int slot, int C, int H, int W, int noise_dim, int tanh_out, const float* blob, size_t n_floats);
int ganrev_forward_G(ganrev_ctx* ctx, const float* noise, int64_t N, float* images);
int ganrev_forward_R(ganrev_ctx* ctx, int slot, const float* images, const uint8_t* mask, int64_t N, float* attrs);
int ganrev_fix_l2(ganrev_ctx* ctx, int slot, const float* images, const uint8_t* mask, int64_t N, float* attrs, float* fixed, double* l2);
int ganrev_l2(ganrev_ctx* ctx, const float* a, const float* b, int64_t N, int px, double* l2);
int ganrev_nearest_l2(ganrev_ctx* ctx, const float* queries, int Q, const float* set, int64_t N, int px, int64_t* ids, double* dist);
int ganrev_anomaly_flags(ganrev_ctx* ctx, const double* l2, int64_t n_calc, int64_t n_show, double quantile, uint8_t* flags, double* thr);
int ganrev_buffer_put(ganrev_ctx* ctx, int which, const void* host, int64_t rows);
int ganrev_buffer_get(ganrev_ctx* ctx, int which, void* host, int64_t row0, int64_t rows);
int ganrev_db_set(ganrev_ctx* ctx, const float* vecs, int64_t N, int d);
int ganrev_cosine(ganrev_ctx* ctx, const float* a, const float* b, int d, float* out);
int ganrev_search_cosine(ganrev_ctx* ctx, const float* queries, int Q, int k, int64_t* ids, float* scores);
int ganrev_search_rows(ganrev_ctx* ctx, const int64_t* rows, int Q, int k, int64_t* ids, float* scores);
int ganrev_kmeans(ganrev_ctx* ctx, int k, int niter, const float* init_centroids, float* centroids, float* total_counts, int32_t* last_labels);
int ganrev_assign_cosine_min(ganrev_ctx* ctx, const float* centroids, int k, int32_t* cluster, float* cosv);
int ganrev_cluster_members(ganrev_ctx* ctx, int k, int m, const float* images, int px, int64_t* member_ids, int32_t* member_counts, float* mean_images);
int ganrev_refine_l2(ganrev_ctx* ctx, int slot, const float* images, const float* z0, int64_t N, int iters, const float* hyper6, float* attrs, float* fixed, double* l2);
int ganrev_train_R_init(ganrev_ctx* ctx, int C, int H, int W, int noise_dim, int tanh_out, int fixer, const float* blob, size_t n_floats);
int ganrev_train_R_step(ganrev_ctx* ctx, const float* noise, int B, const uint8_t* masks, size_t mask_bytes, const float* hyper7, double* loss2);
int ganrev_train_R_state(ganrev_ctx* ctx, int what, float* out, size_t n_floats);
int ganrev_sync(ganrev_ctx* ctx);
int ganrev_set_option(ganrev_ctx* ctx, const char* name, int64_t value);
]]

local lib = ffi.load(os.getenv('GANREV_LIB') or 'ganrev_cuda')   -- libganrev_cuda.so on LD_LIBRARY_PATH
local M = {}

local function check(ctx, rc)
    if rc ~= 0 then error(string.format('ganrev error %d: %s', rc, ffi.string(lib.ganrev_last_error(ctx)))) end
end
local function fptr(t) return t and t:contiguous():data() or nil end   -- FloatTensor:data() -> float*

function M.new(device)
    local out = ffi.new('ganrev_ctx*[1]')
    local rc = lib.ganrev_create(out, device or 0)
    if rc ~= 0 then error('ganrev_create failed (needs an sm_100 GPU; there is no CPU fallback), rc=' .. rc) end
    return ffi.gc(out[0], lib.ganrev_destroy)
end

-- multi-GPU: one Lua state per GPU.  Rank 0 creates the id, the launcher ships the bytes.
function M.unique_id(ctx)
    local buf, len = ffi.new('uint8_t[256]'), ffi.new('size_t[1]')
    check(ctx, lib.ganrev_comm_unique_id(ctx, buf, 256, len))
    return ffi.string(buf, len[0])
end
function M.comm_init(ctx, world, rank, id)
    check(ctx, lib.ganrev_comm_init(ctx, world, rank, id, #id))
end
-- The hand-off as code: one `th apply_r.lua` process per GPU (RANK / WORLD_SIZE in the environment), a path on
-- a file system all of them see.  Rank 0 writes the id to `path .. '.tmp'` and renames it (atomic on POSIX), the
-- others poll for `path`; every rank then joins the communicator.  gan-reverser_b200/dist.py has the same protocol.
function M.comm_init_file(ctx, world, rank, path, timeout_s)
    if world == 1 then return end
    local id
    if rank == 0 then
        id = M.unique_id(ctx)
        local f = assert(io.open(path .. '.tmp', 'wb'))
        f:write(id); f:close()
        assert(os.rename(path .. '.tmp', path))
    else
        local t0 = os.time()
        while true do
            local f = io.open(path, 'rb')
            if f then
                id = f:read('*a'); f:close()
                if #id > 0 then break end
            end
            if os.time() - t0 > (timeout_s or 120) then error('no NCCL unique id at ' .. path) end
            ffi.C.usleep(20000)
        end
    end
    M.comm_init(ctx, world, rank, id)
end

-- Flatten a trained nn.Sequential into the weight blob of include/ganrev.h: every Linear /
-- (cudnn.)SpatialConvolution as weight then bias, every (Spatial)BatchNormalization as
-- gamma, beta, running_mean, running_var -- in module order (models.lua:115-132, 409-451).
function M.flatten(model)
    local parts, n = {}, 0
    local function push(t) t = t:float():contiguous():view(-1); table.insert(parts, t); n = n + t:nElement() end
    for _, m in ipairs(model.modules) do
        local tn = torch.typename(m)
        if tn == 'nn.Linear' or tn:find('SpatialConvolution') then
            push(m.weight); push(m.bias)
        elseif tn:find('BatchNormalization') then
            push(m.weight); push(m.bias); push(m.running_mean)
            -- newer nn keeps running_var, cudnn R3-era nn kept running_std = 1/sqrt(var+eps)
            if m.running_var then push(m.running_var)
            else push(torch.pow(m.running_std:float(), -2):add(-(m.eps or 1e-5))) end
        end
    end
    local blob, o = torch.FloatTensor(n), 1
    for _, t in ipairs(parts) do blob:narrow(1, o, t:nElement()):copy(t); o = o + t:nElement() end
    return blob
end

-- Weight blobs without nn / cudnn -----------------------------------------------------------
-- Layout of include/ganrev.h ("Weight blob"), as {kind, n_out, fan_in} records in models.lua module order.
local function g_layout(C, H, W, nd)
    local F = 512 * (H / 4) * (W / 4)
    return {{'w', F, nd}, {'bn', F}, {'w', 256, 512 * 9}, {'bn', 256}, {'w', 128, 256 * 9}, {'bn', 128}, {'w', C, 128 * 9}}
end
local function r_layout(C, H, W, nd)
    local F = 128 * (H / 4) * (W / 4)
    return {{'w', 64, C * 9}, {'bn', 64}, {'w', 64, 64 * 9}, {'bn', 64}, {'w', 64, 64 * 9}, {'bn', 64}, {'w', 128, 64 * 9}, {'bn', 128},
            {'w', 128, 128 * 9}, {'bn', 128}, {'w', 128, 128 * 9}, {'bn', 128}, {'w', 512, F}, {'bn', 512}, {'w', nd, 512}}
end
-- Random init = what models.lua + w_init(net, 'heuristic') leave behind (weight-init.lua:14-16, 52-73): weights
-- U(+-1/sqrt(fan_in)), every bias (BN beta included) zero, BN gamma U(0,1), running mean 0 / var 1.  Drawn from
-- torch's global generator, so torch.manualSeed(OPT.seed) (apply_r.lua:35) makes it reproducible.
local function init_blob(layout)
    local n = 0
    for _, l in ipairs(layout) do n = n + (l[1] == 'w' and l[2] * l[3] + l[2] or 4 * l[2]) end
    local blob, o = torch.FloatTensor(n):zero(), 1
    for _, l in ipairs(layout) do
        if l[1] == 'w' then
            local bound = 1 / math.sqrt(l[3])
            blob:narrow(1, o, l[2] * l[3]):uniform(-bound, bound); o = o + l[2] * l[3] + l[2]      -- bias stays zero
        else
            blob:narrow(1, o, l[2]):uniform(0, 1)                                                -- gamma
            blob:narrow(1, o + 3 * l[2], l[2]):fill(1); o = o + 4 * l[2]                          -- running_var
        end
    end
    return blob
end
function M.init_blob_G(dimensions, noiseDim) return init_blob(g_layout(dimensions[1], dimensions[2], dimensions[3], noiseDim)) end
function M.init_blob_R(dimensions, noiseDim) return init_blob(r_layout(dimensions[1], dimensions[2], dimensions[3], noiseDim)) end
-- A trained checkpoint converted offline by `python tools/net2blob.py logs/adversarial.net` (Torch7 .net -> raw float32
-- blob + a .json with the geometry): the Lua process then needs neither nn nor cudnn to deserialise it.
function M.read_blob(path)
    return torch.FloatTensor(torch.FloatStorage(path))
end

-- MODELS.create_G(dimensions, noiseDim, cuda)   models.lua:201-203: random-init G3 living in the library
function M.create_G(ctx, dimensions, noiseDim, blob)
    return M.wrap_G(ctx, blob or M.init_blob_G(dimensions, noiseDim), dimensions, noiseDim)
end
-- MODELS.create_R(dimensions, noiseDim, noiseMethod, fixer, cuda)   models.lua:385-387
function M.create_R(ctx, dimensions, noiseDim, noiseMethod, fixer, blob)
    return M.wrap_R(ctx, blob or M.init_blob_R(dimensions, noiseDim), fixer and 1 or 0, dimensions, noiseDim, noiseMethod, fixer)
end

-- Object with the nn.Module protocol apply_r.lua uses (:forward, :evaluate, :training, :float) over a trained
-- nn.Sequential (flattened here) or a ready weight blob (a torch.FloatTensor).
function M.wrap_G(ctx, model, dimensions, noiseDim)
    local blob = torch.isTensor(model) and model:float():contiguous() or M.flatten(model)
    check(ctx, lib.ganrev_load_G(ctx, dimensions[1], dimensions[2], dimensions[3], noiseDim, blob:data(), blob:nElement()))
    local G = {ctx = ctx, dimensions = dimensions, noiseDim = noiseDim}
    function G:forward(noise)                                  -- utils/nn_utils.lua:5-33 batches; the library chunks internally
        noise = noise:float():contiguous()
        if noise:dim() == 1 then noise = noise:view(1, -1) end
        local N = noise:size(1)
        local images = torch.FloatTensor(N, dimensions[1], dimensions[2], dimensions[3])
        check(ctx, lib.ganrev_forward_G(ctx, noise:data(), N, images:data()))
        self.output = images
        return images
    end
    function G:evaluate() return self end
    function G:training() error('libganrev_cuda implements inference only') end
    function G:float() error('no CPU fallback: the apply_r path runs on the B200 only') end
    function G:cuda() return self end
    return G
end

-- MODELS.create_R(dimensions, noiseDim, noiseMethod, fixer, cuda) replacement.  slot 0 = R,
-- slot 1 = R_fixer.  The fixer's always-on input Dropout(0.5) (models.lua:399-406) is drawn
-- here with torch.bernoulli and passed down as an explicit mask (x*mask, no rescale).
function M.wrap_R(ctx, model, slot, dimensions, noiseDim, noiseMethod, fixer)
    assert(noiseMethod == 'normal' or noiseMethod == 'uniform')          -- models.lua:390
    local blob = torch.isTensor(model) and model:float():contiguous() or M.flatten(model)
    check(ctx, lib.ganrev_load_R(ctx, slot, dimensions[1], dimensions[2], dimensions[3], noiseDim,
                                 noiseMethod ~= 'normal' and 1 or 0, blob:data(), blob:nElement()))
    local R = {ctx = ctx, slot = slot, fixer = fixer, noiseDim = noiseDim}
    function R:forward(images, mask)
        images = images:float():contiguous()
        if images:dim() == 3 then images = images:view(1, images:size(1), images:size(2), images:size(3)) end
        local N = images:size(1)
        if self.fixer and mask == nil then
            mask = torch.ByteTensor(images:size()):bernoulli(0.5)
        end
        local attrs = torch.FloatTensor(N, noiseDim)
        check(ctx, lib.ganrev_forward_R(ctx, slot, images:data(), mask and mask:contiguous():data() or nil, N, attrs:data()))
        self.output = attrs
        return attrs
    end
    function R:evaluate() return self end
    function R:training() error('libganrev_cuda implements inference only') end
    function R:float() error('no CPU fallback: the apply_r path runs on the B200 only') end
    function R:cuda() return self end
    return R
end

-- cosineSimilarity(v1, v2)  apply_r.lua:396-400
function M.cosineSimilarity(ctx, v1, v2)
    local out = ffi.new('float[1]')
    v1, v2 = v1:float():contiguous(), v2:float():contiguous()
    check(ctx, lib.ganrev_cosine(ctx, v1:data(), v2:data(), v1:nElement(), out))
    return tonumber(out[0])
end

-- unsup.kmeans(x, k, niter)  apply_r.lua:198 -> centroids, counts.  The N(0,1) row-normalised
-- initial centroids unsup draws internally are drawn here (same torch RNG stream position).
function M.kmeans(ctx, x, k, niter, init)
    x = x:float():contiguous()
    local N, d = x:size(1), x:size(2)
    if not init then
        init = torch.FloatTensor(k, d):normal()
        for i = 1, k do init[i]:div(init[i]:norm()) end
    end
    check(ctx, lib.ganrev_db_set(ctx, x:data(), N, d))
    local cen, counts = torch.FloatTensor(k, d), torch.FloatTensor(k)
    check(ctx, lib.ganrev_kmeans(ctx, k, niter, init:contiguous():data(), cen:data(), counts:data(), nil))
    return cen, counts
end

-- createClusterImages inner loops  apply_r.lua:206-243.  Returns 1-based img2cluster, the
-- per-cluster member lists (1-based, sorted by cosine descending) and the mean faces.
function M.cluster(ctx, attributes, centroids, images, nbMaxPerCluster)
    attributes, images = attributes:float():contiguous(), images:float():contiguous()
    local N, k = attributes:size(1), centroids:size(1)
    check(ctx, lib.ganrev_db_set(ctx, attributes:data(), N, attributes:size(2)))
    local cl, cv = torch.IntTensor(N), torch.FloatTensor(N)
    check(ctx, lib.ganrev_assign_cosine_min(ctx, centroids:float():contiguous():data(), k, cl:data(), cv:data()))
    local px = images:nElement() / N
    local ids, cnt = torch.LongTensor(k, nbMaxPerCluster), torch.IntTensor(k)
    local mean = torch.FloatTensor(k, px)
    check(ctx, lib.ganrev_cluster_members(ctx, k, nbMaxPerCluster, images:data(), px, ids:data(), cnt:data(), mean:data()))
    return cl:add(1), cv, ids:add(1), cnt, mean
end

-- createSimilaritySearchImages inner loops  apply_r.lua:267-282: ids (1-based) and scores of the
-- k most similar database rows for each query row.
function M.search(ctx, db, queries, k)
    db, queries = db:float():contiguous(), queries:float():contiguous()
    check(ctx, lib.ganrev_db_set(ctx, db:data(), db:size(1), db:size(2)))
    local Q = queries:size(1)
    local ids, scores = torch.LongTensor(Q, k), torch.FloatTensor(Q, k)
    check(ctx, lib.ganrev_search_cosine(ctx, queries:data(), Q, k, ids:data(), scores:data()))
    return ids:add(1), scores
end

-- the same with the needles given as (1-based) rows of db itself, apply_r.lua:268
function M.search_rows(ctx, db, needle_rows, k)
    db = db:float():contiguous()
    check(ctx, lib.ganrev_db_set(ctx, db:data(), db:size(1), db:size(2)))
    local Q = needle_rows:size(1)
    local rows0 = needle_rows:long():add(-1):contiguous()
    local ids, scores = torch.LongTensor(Q, k), torch.FloatTensor(Q, k)
    check(ctx, lib.ganrev_search_rows(ctx, rows0:data(), Q, k, ids:data(), scores:data()))
    return ids:add(1), scores
end

-- detectAnomalies  apply_r.lua:355-378: fixed = G(attributesFixer); dist = torch.dist per image;
-- flags = (1 - dist) <= sorted[floor(n*threshold)]
function M.anomalies(ctx, images, fixed, nbImagesCalculations, nbImagesShow, threshold)
    images, fixed = images:float():contiguous(), fixed:float():contiguous()
    local n = nbImagesCalculations
    local px = images:nElement() / images:size(1)
    local l2 = torch.DoubleTensor(n)
    check(ctx, lib.ganrev_l2(ctx, images:data(), fixed:data(), n, px, l2:data()))
    local flags, thr = torch.ByteTensor(nbImagesShow), ffi.new('double[1]')
    check(ctx, lib.ganrev_anomaly_flags(ctx, l2:data(), n, nbImagesShow, threshold, flags:data(), thr))
    return flags, l2:mul(-1):add(1), tonumber(thr[0])
end

-- New work (the reference stops at R's single pass, apply_r.lua:152-153): refine recovered vectors by gradient descent through G.
-- images = N x C x H x W, attributes = N x noiseDim (R's or R_fixer's output, the starting point), nbIterations Adam steps on
-- ||G(z) - x||^2 + prior ||z||^2 per image; opt = {lr, beta1, beta2, eps, prior, zclamp} (defaults 0.01, 0.9, 0.999, 1e-8, 0, 0 = no
-- clamp).  slot = which ATTRS buffer keeps the result (default 1, the fixer's).  Returns refined attributes, G(refined), distances.
function M.refine_l2(ctx, images, attributes, nbIterations, opt, slot)
    opt = opt or {}
    images, attributes = images:float():contiguous(), attributes:float():contiguous()
    local N = images:size(1)
    local hyper = torch.FloatTensor({opt.lr or 0.01, opt.beta1 or 0.9, opt.beta2 or 0.999, opt.eps or 1e-8, opt.prior or 0, opt.zclamp or 0})
    local refined, fixed, l2 = torch.FloatTensor(N, attributes:size(2)), torch.FloatTensor(images:size()), torch.DoubleTensor(N)
    check(ctx, lib.ganrev_refine_l2(ctx, slot or 1, images:data(), attributes:data(), N, nbIterations, hyper:data(),
                                    refined:data(), fixed:data(), l2:data()))
    return refined, fixed, l2
end

-- findClosestNeighboursOf  sample.lua:128-148: images = list of image tensors, trainingSet = N x C x H x W tensor.
-- Returns the same list of {image, closest training image, distance}.
function M.findClosestNeighboursOf(ctx, images, trainingSet)
    local Q = #images
    if Q == 0 then return {} end
    local q = torch.FloatTensor(Q, images[1]:nElement())
    for i = 1, Q do q[i]:copy(images[i]:float():view(-1)) end
    local ts = trainingSet:float():contiguous()
    local N, px = ts:size(1), ts:nElement() / ts:size(1)
    local ids, dist = torch.LongTensor(Q), torch.DoubleTensor(Q)
    check(ctx, lib.ganrev_nearest_l2(ctx, q:data(), Q, ts:data(), N, px, ids:data(), dist:data()))
    local result = {}
    for i = 1, Q do
        table.insert(result, {images[i], ts[ids[i] + 1]:clone(), dist[i]})
    end
    return result
end

-- train_r.lua:129-170.  trainer = ganrev.train_R(ctx, dimensions, noiseDim, noiseMethod, fixer, blob): the optimiser state (Adam's
-- m / v, step count) lives in the context; G must be loaded (train_r.lua:96-98).  trainer.step(noise, masks, hyper) replaces
--   optim.adam(fevalR, PARAMETERS_R, OPTSTATE.adam.R)   train_r.lua:165
-- noise = NN_UTILS.createNoiseInputs(OPT.batchSize); masks = list of ByteTensors in module order (include/ganrev.h), drawn by the
-- caller with torch.bernoulli so Torch's generator keeps owning the randomness; hyper = {learningRate, beta1, beta2, epsilon,
-- R_L1, R_L2, R_clamp} (defaults: optim.adam's + train_r.lua:22-24).  Returns the criterion's loss and feval's f (with penalties).
function M.train_R(ctx, dimensions, noiseDim, noiseMethod, fixer, blob)
    blob = (blob or M.init_blob_R(dimensions, noiseDim)):float():contiguous()
    check(ctx, lib.ganrev_train_R_init(ctx, dimensions[1], dimensions[2], dimensions[3], noiseDim,
                                       noiseMethod ~= 'normal' and 1 or 0, fixer and 1 or 0, blob:data(), blob:nElement()))
    local n_floats = blob:nElement()
    local T = {}
    function T.step(noise, masks, hyper)
        local z = noise:float():contiguous()
        local total = 0
        for _, m in ipairs(masks) do total = total + m:nElement() end
        local mk = torch.ByteTensor(total)
        local at = 1
        for _, m in ipairs(masks) do mk:narrow(1, at, m:nElement()):copy(m:byte():view(-1)); at = at + m:nElement() end
        local hy = torch.FloatTensor(hyper or {1e-3, 0.9, 0.999, 1e-8, 0, 1e-4, 1})
        local out = ffi.new('double[2]')
        check(ctx, lib.ganrev_train_R_step(ctx, z:data(), z:size(1), mk:data(), total, hy:data(), out))
        return tonumber(out[0]), tonumber(out[1])
    end
    -- what: 0 parameters + running statistics (the blob create_R / ganrev_load_R take, what train_r.lua:228-235 saves),
    -- 1 last gradients, 2 / 3 Adam's m / v
    function T.state(what)
        local out = torch.FloatTensor(n_floats)
        check(ctx, lib.ganrev_train_R_state(ctx, what or 0, out:data(), n_floats))
        return out
    end
    return T
end

return M
